#!/usr/bin/env python
"""Generate the golden fixtures of tests/golden/ by running THE REFERENCE'S OWN CUDA KERNELS (oracle/_ref, built from a checkout
of the reference by oracle/build_ref.py for sm_100a) on seeded inputs.  Run on a B200:

    python tests/golden/make_golden.py OUTDIR      # then copy OUTDIR/*.npz to tests/golden/

Inputs are regenerated from seeds by the tests (tests/_golden_inputs.py); only outputs (and tiny inputs) are stored, so the
fixtures stay small.  The reference has no golden vectors or tests of its own (SURVEY.md section 4); these files are what
pins the CPU oracle (tests/test_oracle_cpu.py compares oracle/ntx_oracle.c against them without any GPU).

tests/golden/reference_outputs.npz, what the GPU tests compare with the reference's kernels, is written by those tests themselves
(tests/_util.py: reference_output), on a B200 with oracle/_ref built:

    NTX_RECORD_REFERENCE=$PWD/tests/golden/reference_outputs.npz python -m pytest -m gpu \
        tests/test_gpu_grid.py tests/test_gpu_mlp.py tests/test_gpu_training.py tests/test_gpu_field.py tests/test_gpu_sh.py tests/test_gpu_raymarching.py
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from _golden_inputs import GRID_CASES, MLP_CASES, grid_case_inputs, mlp_case_inputs, scene_inputs, sh_inputs  # noqa: E402
from _util import _digest, ref  # noqa: E402

DEV = "cuda"
SAMPLE = 512


def shrink_grid(out, name):
    """keep grid.npz small: the outputs as a digest of the whole array plus a fixed seeded sample of its elements, the table and
    input gradients as a seeded sample of rows plus the largest magnitude of the whole"""
    rng = np.random.default_rng(0)
    for k in ("_out_LBC", "_dy_dx"):
        a = out.pop(name + k).reshape(-1)
        a = a.view({2: np.uint16, 4: np.uint32}[a.itemsize])          # compared bit for bit
        idx = np.sort(rng.choice(a.size, SAMPLE, replace=False))
        out[name + k + ":rows"], out[name + k + ":sample"], out[name + k + ":digest"] = idx.astype(np.int32), a[idx], _digest(a)
    rows, vals = out.pop(name + "_grad_rows"), out.pop(name + "_grad_vals")
    sel = np.sort(rng.choice(len(rows), min(SAMPLE, len(rows)), replace=False))
    out[name + "_grad_rows"], out[name + "_grad_vals"] = rows[sel].astype(np.int32), vals[sel]
    out[name + "_grad_vals_absmax"] = np.abs(vals.astype(np.float64)).max()
    gi = out.pop(name + "_grad_inputs")
    sel = np.sort(rng.choice(len(gi), min(SAMPLE, len(gi)), replace=False))
    out[name + "_grad_inputs:rows"], out[name + "_grad_inputs:sample"] = sel.astype(np.int32), gi[sel]
    out[name + "_grad_inputs_absmax"] = np.abs(gi.astype(np.float64)).max()


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def main(outdir):
    os.makedirs(outdir, exist_ok=True)
    g, f, s, r = ref("gridencoder"), ref("ffmlp"), ref("shencoder"), ref("raymarching")

    # ---- the device's per-level scales (exp2f is an approximate instruction on the GPU) ---------------------------
    import nerf_texture_b200
    from nerf_texture_b200 import _lib as L
    out = {}
    for name, case in GRID_CASES.items():
        x, emb, offsets, pls, cfg = grid_case_inputs(case)
        nlev = offsets.shape[0] - 1
        sc = torch.empty(nlev, device=DEV)
        L.call("ntx_grid_level_scales", float(np.log2(pls)), cfg["base_resolution"], nlev, sc.data_ptr(), L.stream())
        B, D = x.shape
        C = emb.shape[1]
        xt, et, ot = T(x), T(emb), T(offsets)
        o = torch.empty(nlev, B, C, dtype=et.dtype, device=DEV)
        dy = torch.empty(B, nlev * D * C, dtype=et.dtype, device=DEV)
        g.grid_encode_forward(xt, et, ot, o, B, D, C, nlev, float(np.log2(pls)), cfg["base_resolution"], True, dy, case["gridtype"], cfg["align_corners"])
        grad = T(np.random.default_rng(case["seed"] + 100).standard_normal((nlev, B, C)).astype(emb.dtype))
        ge = torch.zeros_like(et)
        gi = torch.zeros(B, D, dtype=et.dtype, device=DEV)
        g.grid_encode_backward(grad, xt, et, ot, ge, B, D, C, nlev, float(np.log2(pls)), cfg["base_resolution"], True, dy, gi, case["gridtype"], cfg["align_corners"])
        torch.cuda.synchronize()
        out[name + "_scales"] = sc.cpu().numpy()
        out[name + "_out_LBC"] = o.cpu().numpy()
        out[name + "_dy_dx"] = dy.cpu().numpy()
        nz = torch.nonzero(ge.float().abs().sum(1)).flatten().cpu().numpy()[:4096]      # sparse sample of the table gradient
        out[name + "_grad_rows"] = nz.astype(np.int64)
        out[name + "_grad_vals"] = ge[torch.from_numpy(nz).to(DEV)].cpu().numpy()
        out[name + "_grad_inputs"] = gi.cpu().numpy()
        shrink_grid(out, name)
    np.savez_compressed(os.path.join(outdir, "grid.npz"), **out)

    out = {}
    for name, case in MLP_CASES.items():
        x, w = mlp_case_inputs(case)
        B = x.shape[0]
        f.allocate_splitk(case["layers"] + 1)
        o = torch.empty(B, 16, dtype=torch.half, device=DEV)
        buf = torch.empty(B, case["hidden"], dtype=torch.half, device=DEV)
        f.ffmlp_inference(T(x), T(w), B, case["in_dim"], 16, case["hidden"], case["layers"], 0, 6, buf, o)
        fb = torch.empty(case["layers"], B, case["hidden"], dtype=torch.half, device=DEV)
        o2 = torch.empty(B, 16, dtype=torch.half, device=DEV)
        f.ffmlp_forward(T(x), T(w), B, case["in_dim"], 16, case["hidden"], case["layers"], 0, 6, fb, o2)
        torch.cuda.synchronize()
        out[name + "_out"] = o.cpu().numpy()
        out[name + "_fwd_last"] = fb[-1].cpu().numpy()
    np.savez_compressed(os.path.join(outdir, "ffmlp.npz"), **out)

    out = {}
    for deg in (1, 2, 4, 6, 8):
        d = sh_inputs(deg)
        B = d.shape[0]
        o = torch.empty(B, deg * deg, device=DEV)
        dy = torch.empty(B, 3 * deg * deg, device=DEV)
        s.sh_encode_forward(T(d), o, B, 3, deg, True, dy)
        torch.cuda.synchronize()
        out["deg%d_out" % deg] = o.cpu().numpy()
        out["deg%d_dy_dx" % deg] = dy.cpu().numpy()
    np.savez_compressed(os.path.join(outdir, "sh.npz"), **out)

    out = {}
    for name in ("c1", "c2"):
        sc = scene_inputs(name)
        o, d, bits, aabb = T(sc["rays_o"]), T(sc["rays_d"]), T(sc["bits"]), T(sc["aabb"])
        N = sc["rays_o"].shape[0]
        nears, fars = torch.empty(N, device=DEV), torch.empty(N, device=DEV)
        r.near_far_from_aabb(o, d, aabb, N, 0.2, nears, fars)
        M = N * sc["max_steps"]
        xyzs, dirs, deltas = torch.zeros(M, 3, device=DEV), torch.zeros(M, 3, device=DEV), torch.zeros(M, 2, device=DEV)
        rays = torch.empty(N, 3, dtype=torch.int32, device=DEV)
        cnt = torch.zeros(2, dtype=torch.int32, device=DEV)
        r.march_rays_train(o, d, bits, sc["bound"], sc["dt_gamma"], sc["max_steps"], N, sc["cascade"], sc["H"], M, nears, fars, xyzs, dirs, deltas, rays, cnt, sc["perturb"])
        torch.cuda.synchronize()
        rays_np = rays.cpu().numpy()
        order = np.argsort(rays_np[:, 0], kind="stable")     # the reference's row order is arbitrary (atomics): store sorted by ray id
        m = int(cnt[0].item())
        rng = np.random.default_rng(7)
        sig = (rng.random(m + 128).astype(np.float32) * 20)
        rgb = rng.random((m + 128, 3)).astype(np.float32)
        ws, dp, im = torch.empty(N, device=DEV), torch.empty(N, device=DEV), torch.empty(N, 3, device=DEV)
        r.composite_rays_train_forward(T(sig), T(rgb), deltas[:m + 128].contiguous(), rays, m + 128, N, ws, dp, im)
        torch.cuda.synchronize()
        out[name + "_nears"], out[name + "_fars"] = nears.cpu().numpy(), fars.cpu().numpy()
        out[name + "_counter"] = cnt.cpu().numpy()
        out[name + "_ray_counts"] = rays_np[order][:, 2]
        # per-ray samples in ray order (what an ordered allocation produces)
        xs, ds = xyzs.cpu().numpy(), deltas.cpu().numpy()
        segs_x = [xs[a:a + c] for a, c in zip(rays_np[order][:, 1], rays_np[order][:, 2])]
        segs_d = [ds[a:a + c] for a, c in zip(rays_np[order][:, 1], rays_np[order][:, 2])]
        out[name + "_xyzs_ordered"] = np.concatenate(segs_x) if m else np.zeros((0, 3), np.float32)
        out[name + "_deltas_ordered"] = np.concatenate(segs_d) if m else np.zeros((0, 2), np.float32)
        out[name + "_ws"], out[name + "_depth"], out[name + "_image"] = ws.cpu().numpy(), dp.cpu().numpy(), im.cpu().numpy()
        out[name + "_comp_ray_order"] = rays_np[:, 0]         # which image row each reference ray row wrote (needed to re-index sig/rgb)
        out[name + "_comp_offsets"] = rays_np[:, 1]
        # one inference-loop iteration: march_rays (n_step 4) + composite_rays + compact_rays
        alive = torch.arange(N, dtype=torch.int32, device=DEV)
        tt = nears.clone()
        n_step = 4
        Mi = N * n_step + 128 - (N * n_step) % 128
        ix, idr, idl = torch.zeros(Mi, 3, device=DEV), torch.zeros(Mi, 3, device=DEV), torch.zeros(Mi, 2, device=DEV)
        r.march_rays(N, n_step, alive, tt, o, d, sc["bound"], sc["dt_gamma"], sc["max_steps"], sc["cascade"], sc["H"], bits, nears, fars, ix, idr, idl, sc["perturb"])
        sig2 = T(rng.random(Mi).astype(np.float32) * 200)
        rgb2 = T(rng.random((Mi, 3)).astype(np.float32))
        ws2, dp2, im2 = torch.zeros(N, device=DEV), torch.zeros(N, device=DEV), torch.zeros(N, 3, device=DEV)
        r.composite_rays(N, n_step, alive, tt, sig2, rgb2, idl, ws2, dp2, im2)
        alive2, t2 = torch.zeros_like(alive), torch.zeros_like(tt)
        c2 = torch.zeros(1, dtype=torch.int32, device=DEV)
        r.compact_rays(N, alive2, alive, t2, tt, c2)
        torch.cuda.synchronize()
        k = int(c2.item())
        a2, t2n = alive2[:k].cpu().numpy(), t2[:k].cpu().numpy()
        o2 = np.argsort(a2, kind="stable")
        out[name + "_inf_xyzs"], out[name + "_inf_deltas"] = ix.cpu().numpy(), idl.cpu().numpy()
        out[name + "_inf_t_after"] = tt.cpu().numpy()
        out[name + "_inf_ws"], out[name + "_inf_image"], out[name + "_inf_depth"] = ws2.cpu().numpy(), im2.cpu().numpy(), dp2.cpu().numpy()
        out[name + "_inf_alive_sorted"], out[name + "_inf_t_sorted"] = a2[o2], t2n[o2]
    np.savez_compressed(os.path.join(outdir, "raymarching.npz"), **out)
    for fn in sorted(os.listdir(outdir)):
        print(fn, os.path.getsize(os.path.join(outdir, fn)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE))
