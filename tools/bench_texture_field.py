#!/usr/bin/env python
"""Fused texture-field density (ntx_texture_field_density) against the same computation composed from the in-tree drop-ins:

    python tools/bench_texture_field.py [--lat 340] [--iters 10]

Two workloads on the 230 K-triangle bumpy sphere of tools/bench_mesh.py, bound 1, cfgT texture grid, the tinycudann shim's sigma_net
(41 -> 32 -> 16), h_threshold 0.1, under fp16 autocast without gradients (how update_extra_state calls NeRFNetwork.density):
  (a) `shell`: 2^20 samples of 8192 camera-like rays x 128 steps through 0.45 <= |x| <= 0.95, in ray order (bench_mesh.py's generator);
  (b) `grid`: the 128^3 cell centres of a full density-grid update of cascade 0 (renderer.py:585-600: 2 * coords / (H - 1) - 1, scaled
      by bound - half_grid_size), in one call — the renderer's chunk S = 128 covers the whole 128^3 grid.
Arms: `composed` = Mesh.project -> GridEncoder -> frequency encoding -> tinycudann.Network -> exp / where; `fused` = texture.density.
Both visit batches of mesh.SORT_MIN samples or more in Morton order.  CUDA events, 3 warm-up calls, a 256 MB write between timed calls
flushes L2, the two arms alternate, median of --iters.  The outputs of both arms are compared bit for bit at the timed size.  Prints
`RESULT {json}` with the GPU's name and power limit.  Reads nothing outside this repository."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _gpu():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in q.stdout.strip().split(",")]
        return name, power
    except Exception as e:                                    # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(e).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lat", type=int, default=340)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--log2-samples", type=int, default=20)
    args = ap.parse_args()
    import numpy as np
    import torch
    import _util as U
    import nerf_texture_b200
    nerf_texture_b200.install()
    from nerf_texture_b200 import texture
    from test_gpu_texture_field import Field, Model, Projector
    assert torch.cuda.is_available(), "this benchmark needs a GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)

    v, f, vn = U.bumpy_sphere(args.lat, args.lat)
    model = Model(Field(Projector(v, f, vn)))

    # (a) shell samples in ray order (tools/bench_mesh.py)
    N = 1 << args.log2_samples
    steps = 128
    rays = N // steps
    g = torch.Generator(device="cpu").manual_seed(0)
    o = torch.nn.functional.normalize(torch.randn(rays, 3, generator=g), dim=-1) * 1.5
    tgt = torch.nn.functional.normalize(torch.randn(rays, 3, generator=g), dim=-1) * 0.6
    d = torch.nn.functional.normalize(tgt - o, dim=-1)
    ts = torch.linspace(0.4, 2.4, steps)
    x = (o[:, None] + ts[None, :, None] * d[:, None]).reshape(-1, 3)
    rad = x.norm(dim=-1)
    shell = torch.where(((rad < 0.45) | (rad > 0.95))[:, None], x / rad[:, None] * rad.clamp(0.45, 0.95)[:, None], x).contiguous().to(dev)
    # (b) cell centres of cascade 0 of a 128^3 density grid, bound 1 (renderer.py:585-598, no jitter)
    H, bound = 128, 1.0
    c = torch.arange(H, dtype=torch.int32, device=dev)
    X, Y, Z = torch.meshgrid(c, c, c, indexing="ij")
    coords = torch.stack([X.reshape(-1), Y.reshape(-1), Z.reshape(-1)], -1)
    hgs = bound / H
    cells = ((2 * coords.float() / (H - 1) - 1) * (bound - hgs)).contiguous()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    arms = {"composed": lambda q: model.density(q), "fused": lambda q: texture.density(model, q)}
    result = {}
    name, power = _gpu()
    with torch.no_grad(), torch.autocast("cuda", torch.float16):
        for wl, q in (("shell", shell), ("grid", cells)):
            outs = {}
            for arm, fn in arms.items():
                for _ in range(3):
                    outs[arm] = fn(q)
            torch.cuda.synchronize()
            assert model.calls > 0
            same = (torch.equal(outs["fused"]["sigma"].view(torch.int32), outs["composed"]["sigma"].view(torch.int32))
                    and torch.equal(outs["fused"]["geo_feat"].view(torch.int16), outs["composed"]["geo_feat"].view(torch.int16)))
            ms = {a: [] for a in arms}
            for _ in range(args.iters):
                for arm, fn in arms.items():
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn(q)
                    e1.record()
                    torch.cuda.synchronize()
                    ms[arm].append(e0.elapsed_time(e1))
            med = {a: float(np.median(t)) for a, t in ms.items()}
            result[wl] = {"samples": int(q.shape[0]), "composed_ms": med["composed"], "fused_ms": med["fused"],
                          "fused_over_composed": med["fused"] / med["composed"], "outputs_equal": bool(same),
                          "in_shell": float((outs["fused"]["sigma"] > 0).float().mean().item()),
                          "composed_ms_all": [round(t, 4) for t in ms["composed"]], "fused_ms_all": [round(t, 4) for t in ms["fused"]]}
            print("%-6s N=%-8d composed %.3f ms  fused %.3f ms  fused/composed %.3f  outputs equal: %s" % (
                wl, q.shape[0], med["composed"], med["fused"], med["fused"] / med["composed"], same), flush=True)
    result.update({"gpu": name, "power_limit": power, "mesh_triangles": int(len(f)), "iters": args.iters})
    print("RESULT " + json.dumps(result))


if __name__ == "__main__":
    main()
