#!/usr/bin/env python
"""bench.py — ray-samples/sec of the per-ray-sample hot path (march -> hash-grid -> fused MLPs -> composite) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one 1024x1024 frame of BASELINE config 3 (random-weight network_ff field, ball occupancy, bound 1, dt_gamma 0,
max_steps 1024) rendered through the libntx C ABI; with N > 1 the frame's rays are sharded over the ranks in interleaved
tiles and the result is all-gathered (config 4, strong scaling).  `value` = non-sentinel samples of the frame / device
time (CUDA events, max over ranks, inputs resident in HBM); `e2e` = the same with rays coming from pinned host memory and
the image read back every step.  `roofline` is for the dominant kernel (the fused field kernel: hash-grid gather + both
MLPs), measured live with CUDA events around every launch of one extra frame.  `cfg2` reports BASELINE config 2 (2^20
random and ray-coherent samples through the fused field kernel and through the stand-alone grid encoder).
`cpu_baseline` / `--impl reference`: the reference has no CPU implementation of this path (SURVEY F1), so the CPU arm is
the oracle port (oracle/ntx_oracle.c, OpenMP over all host cores) rendering a strided sub-sample of the same frame.
`--dump-outputs DIR` writes the frame the last timed step returned (image, depth, weights_sum) as DIR/<name>.npy in float32; the
scene is seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ray-samples/sec (encoder+MLP+composite)"
UNIT = "samples/s"
IMG = 1024
FIELD_BYTES_PER_SAMPLE = 12 + 12 + 4 + 512 + 4 + 12   # xyz, dir, delta | 16 levels x 8 corners x 2 x fp16 | sigma, rgb  (DESIGN.md)
GRID_BYTES_PER_SAMPLE = 12 + 512 + 64                 # SURVEY.md 8d: stand-alone encoder, fp16 table


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """samples nvidia-smi SM clocks + throttle reasons while the timed region runs"""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        # NVML from a thread (a sample every ~5 ms: a timed region of ten 8 ms frames gets ~16 of them); nvidia-smi -lms as fallback
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.samples, self.mask, self.running = [], 0, True
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))

            def loop():
                while self.running:
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)))
                        self.mask |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if getattr(self, "nvml", None) is not None:
            self.running = False
            self.thread.join(timeout=1)
            bits = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}
            return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(n for n, b in bits.items() if self.mask & b), "samples": len(self.samples), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_scene(device, seed=0):
    from nerf_texture_b200 import render, scene
    field = render.NGPField.random(device, seed=seed)
    rays_o, rays_d = scene.pinhole_rays(IMG, IMG, device)
    bits = scene.ball_bitfield(1, 128, 1.0, device)
    return field, rays_o, rays_d, bits


def cpu_render_sample(stride=5, steps=1, warmup=0):
    """oracle (CPU) render of every `stride`-th pixel row/column of the same frame; returns samples/s and a description"""
    import numpy as np
    from oracle import oracle as O
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _util import ball_density_grid, pinhole_rays
    o, d = pinhole_rays(IMG, IMG)
    sel = np.zeros((IMG, IMG), bool)
    sel[::stride, ::stride] = True
    o, d = np.ascontiguousarray(o[sel.ravel()]), np.ascontiguousarray(d[sel.ravel()])
    bits = O.packbits(ball_density_grid(1, 128, 1.0), 0.5)
    offs, pls = O.grid_offsets(3, 16, 2, base_resolution=16, log2_hashmap_size=19, desired_resolution=2048, align_corners=True)
    rng = np.random.default_rng(1)
    emb = (rng.random((int(offs[-1]), 2), dtype=np.float32) * 2 - 1).astype(np.float16)
    ws = ((rng.random(64 * (32 + 64 + 16), dtype=np.float32) * 2 - 1) * np.sqrt(3 / 64)).astype(np.float16)
    wc = ((rng.random(64 * (32 + 128 + 16), dtype=np.float32) * 2 - 1) * np.sqrt(3 / 64)).astype(np.float16)
    times, ns = [], 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        _, _, _, ns, _ = O.render_rays(o, d, bits, 1, 128, 1.0, emb, offs, pls, 16, ws, wc)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return ns / dt, dt, ns, O.num_threads(), "oracle port (oracle/ntx_oracle.c, OpenMP): every %dth row/column of the 1024x1024 frame = %d rays, %d samples per step" % (stride, o.shape[0], ns)


def reference_arm(args):
    """`--impl reference`: the CPU port of the reference path on the host cores (the reference itself is CUDA-only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # One OpenMP thread per PHYSICAL core, set before libgomp loads: with the default (one per hardware thread, 128 on the GPU
    # box) the oracle's many short parallel regions ran 10x slower than with 64 threads (measured: 34 K vs 321 K samples/s).
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:
        phys = max(1, (os.cpu_count() or 2) // 2)
    os.environ["OMP_NUM_THREADS"] = str(phys)     # torchrun exports OMP_NUM_THREADS=1 for its workers: override it here
    os.environ.setdefault("OMP_PROC_BIND", "false")
    value, dt, ns, cores, sample = cpu_render_sample(stride=5, steps=max(1, args.steps), warmup=min(1, args.warmup))   # same sub-sample as cpu_baseline
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": "render_1024x1024_network_ff_random_weights (BASELINE config 3), CPU sub-sample", "l2": "n/a (CPU)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ntx", choices=["ntx", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the cfg2 / roofline side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed step returned as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    from nerf_texture_b200 import _lib as L
    from nerf_texture_b200 import render

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    W, K = max(args.warmup, 3), args.steps
    # host side of the rank on the GPU's own NUMA node (pinned staging buffers, frame mailbox, launches); undone for the CPU baseline
    prev_affinity = L.bind_host_thread_to_gpu(local_rank)
    L.lib()
    assert L.lib().ntx_device_ok() == 1, "libntx needs a CC 10.x device"

    field, rays_o, rays_d, bits = build_scene(device)
    N = rays_o.shape[0]
    if world > 1:
        idx = render.shard_indices(N, world, rank).to(device)
        my_o, my_d = rays_o[idx].contiguous(), rays_d[idx].contiguous()
    else:
        my_o, my_d = rays_o, rays_d

    n_max = render._shard_plan(N, world, 1024, device)[1] if world > 1 else None
    # config 4's exchange step: NVLink peer reads fused into the assembly kernel when symmetric memory is available (NTX_EXCHANGE=nccl
    # forces the all-gather), else ONE NCCL all_gather + the assembly kernel
    exchange = render.PeerFrameExchange.create(N, device=device) if (world > 1 and os.environ.get("NTX_EXCHANGE", "peer") != "nccl") else None
    if world > 1:
        flag = torch.tensor([1 if exchange is not None else 0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)                     # all ranks or none
        if int(flag.item()) == 0:
            exchange = None

    def finish(out):
        if world == 1:
            return out
        if exchange is not None:
            res = exchange.assemble(1.0)
            res["iterations"] = out["iterations"]
            return res
        return render.gather_frame(out, N)

    last = {}

    def step_device():
        # this rank's (resident) shard of the frame, rendered straight into its planar send block, + the exchange and the assembly
        # kernel (config 4); one GPU: the frame
        out = render.render_rays(field, my_o, my_d, bits, 1, 128, block_rows=n_max, cache_mip=True, block_out=exchange.block() if exchange is not None else None)
        last["out"] = finish(out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # samples per frame (untimed, counted once: the scene is deterministic)
    cnt = render.render_rays(field, my_o, my_d, bits, 1, 128, count_samples=True)
    n_local = torch.tensor([cnt["n_samples"]], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(n_local)
    samples_per_frame = int(n_local.item())
    iterations = cnt["iterations"]

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)   # > 126 MB L2

    def timed(fn, steps):
        evs = []
        barrier()
        for _ in range(steps):
            flush.zero_()                      # L2 flush between timed iterations (untimed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            evs.append((e0, e1))
        barrier()
        t = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps         # ms per step, max over ranks

    for _ in range(W):
        step_device()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = L.launches
    ms = timed(step_device, K)
    launches = (L.launches - l0) // K
    clocks = sampler.stop() if rank == 0 else None
    value = samples_per_frame / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in last["out"].items():
            if torch.is_tensor(t):
                np.save(os.path.join(args.dump_outputs, name + ".npy"), t.float().cpu().numpy())
    last.clear()

    # ---- end to end: rays from pinned host memory each step, image + depth read back each step --------------------
    h_o, h_d = my_o.cpu().pin_memory(), my_d.cpu().pin_memory()
    d_o, d_d = torch.empty_like(my_o), torch.empty_like(my_d)
    h_img = torch.empty(N, 3, dtype=torch.float32).pin_memory()
    h_dep = torch.empty(N, dtype=torch.float32).pin_memory()

    def step_e2e():
        d_o.copy_(h_o, non_blocking=True); d_d.copy_(h_d, non_blocking=True)
        out = render.render_rays(field, d_o, d_d, bits, 1, 128, block_rows=n_max, cache_mip=True,       # each rank uploads and renders its own shard
                                 block_out=exchange.block() if exchange is not None else None)
        out = finish(out)
        if rank == 0:
            h_img.copy_(out["image"], non_blocking=True); h_dep.copy_(out["depth"], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    step_e2e()
    ms_e2e = timed(step_e2e, max(3, K // 2))
    e2e = {"value": samples_per_frame / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": int(h_o.numel() * 4 * 2 * world), "d2h_bytes_per_step": int(N * 16)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": "render_1024x1024_network_ff_random_weights (BASELINE config 3%s)" % (("; rays sharded in interleaved 1024-ray tiles + " + ("NVLink peer reads fused into the assembly kernel (symmetric memory)" if exchange is not None else "one NCCL all_gather") + ", config 4") if world > 1 else ""),
                   "field": "hashgrid L=16 T=2^19 F=2 fp16 -> FFMLP(32,16,64,2) -> SH4 -> FFMLP(32,3,64,3)", "rays": N, "samples_per_frame": samples_per_frame,
                   "loop_iterations": iterations, "sample_schedule": "n_step = clamp(32N // n_alive, 1, 256) rounded to 4, walk budget %d, rays that cannot reach an occupied cell dropped before the first march (same image as the reference's clamp(N // n_alive, 1, 8): 43 iterations)" % render.WALK_BUDGET,
                   "max_steps": 1024, "dt_gamma": 0, "occupancy": "ball r=0.5, H=128, 1 cascade (its occupancy mip is built once and cached per bit-field version, like the drop-in march_rays)",
                   "l2": "flushed between timed steps (256 MiB memset)", "parallelism": "ray-sharded x%d" % world,
                   "host": "rank thread bound to the GPU's NUMA node (NVML ideal affinity)" if prev_affinity else "no NUMA binding (NVML unavailable)"},
        "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
    }

    # ---- where a rank's time goes at this N (SCALE runs): march / field kernel sums of one frame (CUDA events inside
    #      ntx_render_rays), the rank's whole shard, and the all-gather + assembly — every rank reports, rank 0 prints
    if world > 1:
        flush.zero_()
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        o = render.render_rays(field, my_o, my_d, bits, 1, 128, time_kernels=True, block_rows=n_max, block_out=exchange.block() if exchange is not None else None)
        ev[1].record()
        finish(o)
        ev[2].record()
        torch.cuda.synchronize()
        mine = torch.tensor([o["march_ms"], o["field_ms"], ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), float(o["iterations"])], dtype=torch.float32, device=device)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        line["per_rank_ms"] = [{"rank": r, "march_ms": round(float(v[0]), 3), "field_ms": round(float(v[1]), 3), "shard_ms": round(float(v[2]), 3),
                                "gather_ms": round(float(v[3]), 3), "iterations": int(v[4])} for r, v in enumerate(allr)]

    if rank == 0 and not args.no_extras:
        peaks, peak_src = measured_peaks()
        # ---- roofline of the dominant kernel: every field launch of one frame bracketed by CUDA events -----------------
        # (ntx_render_rays brackets its own march / field launches with CUDA events on the launching stream when asked to:
        #  same code path, schedule and data as the timed step)
        tk = None
        for _ in range(3):
            flush.zero_()
            o = render.render_rays(field, my_o, my_d, bits, 1, 128, count_samples=True, time_kernels=True)
            if tk is None or o["field_ms"] < tk["field_ms"]:
                tk = o
        kt = tk["field_ms"] * 1e-3
        live = tk["n_samples"]
        nlaunch = tk["iterations"]
        achieved = live * FIELD_BYTES_PER_SAMPLE / kt / 1e9
        # DRAM bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum of ALL field-kernel launches of one frame of this build
        # (one ncu pass, tools/gpu/r2_final.sh -> profiles/r02_field_kernel_traffic.json), divided by the launches that did work
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_field_kernel_traffic.json")))
            traffic = int(tj["dram_bytes_all_field_launches_of_one_frame"] / max(nlaunch, 1))
        except Exception:
            pass
        line["roofline"] = {"bound": "hbm", "kernel": "ngp_field_kernel (hash-grid gather + sigma MLP + SH + colour MLP)", "achieved": achieved,
                            "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_src,
                            "algorithmic_bytes_per_launch": live * FIELD_BYTES_PER_SAMPLE / max(nlaunch, 1),
                            "algorithmic_bytes_per_sample": FIELD_BYTES_PER_SAMPLE, "launches": nlaunch, "avg_launch_us": kt / max(nlaunch, 1) * 1e6,
                            "live_samples": live, "kernel_share_of_step": kt * 1e3 / ms, "march_kernel_ms": tk["march_ms"],
                            "msamples_per_s_in_kernel": live / kt / 1e6,
                            "tensor_note": "36864 FLOP/sample on tcgen05: %.1f TFLOP/s achieved inside the kernel" % (live * 36864 / kt / 1e12)}
        # ---- BASELINE config 1: grid_encode forward L=4 T=2^14 F=2 on 4096 random points — the reference has no CPU path (SURVEY F1), so
        #      the "CPU" number is the oracle port on the host cores; the GPU kernel on the same input next to it
        if prev_affinity:
            os.sched_setaffinity(0, prev_affinity)              # CPU legs (cfg1 here, cpu_baseline below) use every host core; the GPU
        line["cfg1"] = bench_cfg1(torch, L, device)             # side measurements that follow are device-timed
        # ---- BASELINE config 2: 2^20 samples through the fused field kernel and the stand-alone encoder ------------
        line["cfg2"] = bench_cfg2(torch, L, field, device, peaks)
        # ---- the reference's own CUDA kernels (rebuilt for sm_100a, oracle/_ref) on the same frame, when the build is present:
        #      context for the headline only — the contract's reference arm (--impl reference) is the CPU oracle
        if world == 1 and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "_ref_raymarching.so")):
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import compare_ref
                line["reference_cuda"] = compare_ref.main(only_frame=True)
            except Exception as e:      # never let the side measurement break the bench line
                line["reference_cuda"] = {"unavailable": repr(e)[:200]}
        # ---- the drop-in path: the reference's UNMODIFIED nerf/renderer.py + nerf/network_ff.py (baseline/_ref/callers) rendering the
        #      same frame through nerf_texture_b200/compat, next to the same files on the reference's own wrappers + CUDA (oracle/_ref)
        if world == 1:
            line["compat"] = run_tool("run_reference_files.py", [["--backend", "ntx", "--size", str(IMG), "--time", "5"],
                                                                 ["--backend", "ref", "--size", str(IMG), "--time", "5"]], ("ntx", "reference_cuda"), "frame_ms")
            # ---- BASELINE config 5: training step (grid + sigma-MLP forward/backward on 2^18 samples) through the operator API
            line["cfg5"] = run_tool("bench_cfg5.py", [["--backend", "ntx"], ["--backend", "ref"]], ("ntx", "reference_cuda"), "step_ms")
            # ---- SURVEY 8 f3, the mesh front end of the texture field: MeshProjector.project on 2^20 samples — one fused kernel vs the
            #      reference's unmodified torch chain on the drop-in frnn / RayTracer packages vs the CPU restatement
            line["mesh"] = run_tool("bench_mesh.py", [[]], ("ntx",), "project_fused_ms").get("ntx")
        if not args.no_cpu_baseline and world == 1:
            if prev_affinity:
                os.sched_setaffinity(0, prev_affinity)          # the CPU arm uses every host core again
            v, dt, ns, cores, sample = cpu_render_sample(stride=5)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "seconds": dt}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_tool(tool, arg_sets, names, key):
    """run tools/<tool> once per argument set in a subprocess (the two operator stacks cannot share a process: both provide
    `gridencoder`, `ffmlp`, ...), collect its RESULT line; speedup = reference / ntx on `key`"""
    out = {}
    for name, extra in zip(names, arg_sets):
        try:
            r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool)] + extra, capture_output=True, text=True, timeout=900)
            res = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
            out[name] = json.loads(res[0][7:]) if res else {"unavailable": (r.stderr or r.stdout)[-300:]}
        except Exception as e:
            out[name] = {"unavailable": repr(e)[:200]}
    if len(names) < 2:
        return out
    a, b = out.get(names[0], {}), out.get(names[1], {})
    if key in a and key in b and a[key] > 0:
        out["speedup_vs_reference_cuda"] = b[key] / a[key]
    return out


def bench_cfg1(torch, L, device):
    import numpy as np
    from oracle import oracle as O
    offs, pls = O.grid_offsets(3, 4, 2, per_level_scale=2, base_resolution=16, log2_hashmap_size=14, align_corners=False)
    rng = np.random.default_rng(1)
    emb = (rng.random((int(offs[-1]), 2), dtype=np.float32) * 2 - 1).astype(np.float32)
    x = np.random.default_rng(0).random((4096, 3), dtype=np.float32)
    ts = []
    for it in range(55):
        t0 = time.perf_counter()
        O.grid_encode(x, emb, offs, pls, 16, gridtype=0, align_corners=False)
        if it >= 5:
            ts.append(time.perf_counter() - t0)
    cpu_us = statistics.median(ts) * 1e6
    xt, et, ot = torch.from_numpy(x).to(device), torch.from_numpy(emb).to(device), torch.from_numpy(np.asarray(offs, np.int32)).to(device)
    out = torch.empty(4096, 8, device=device)
    fn = lambda: L.call("ntx_grid_encode_forward", L.ptr(xt), L.ptr(et), L.ptr(ot), L.ptr(out), 4096, 3, 2, 4, 1.0, 16, 0, None, 0, 0, L.F32, L.LAYOUT_BLC, L.stream())
    for _ in range(5):
        fn()
    evs = []
    for _ in range(50):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    gpu_us = statistics.median(a.elapsed_time(b) for a, b in evs) * 1e3
    return {"cpu_oracle_port_us": cpu_us, "cpu_threads": O.num_threads(), "ntx_gpu_us": gpu_us, "points": 4096,
            "note": "grid_encode forward, L=4 T=2^14 F=2 fp32 table, median of 50; the CPU arm is the oracle port (no reference CPU path exists)"}


def bench_cfg2(torch, L, field, device, peaks):
    import math
    B = 1 << 20
    g = torch.Generator(device="cpu").manual_seed(0)
    x_rand = (torch.rand(B, 3, generator=g) * 2 - 1).to(device)
    d = torch.randn(B, 3, generator=g)
    d = (d / d.norm(dim=1, keepdim=True)).to(device)
    # ray-coherent variant: 4096 rays x 256 steps of dt_min through the unit cube
    o = (torch.rand(4096, 1, 3, generator=g) * 0.6 - 0.3)
    dd = torch.randn(4096, 1, 3, generator=g); dd = dd / dd.norm(dim=-1, keepdim=True)
    t = (torch.arange(256).float() * (2 * math.sqrt(3) / 1024)).view(1, 256, 1)
    x_coh = (o + dd * t).clamp(-1, 1).reshape(-1, 3).contiguous().to(device)
    d_coh = dd.expand(4096, 256, 3).reshape(-1, 3).contiguous().to(device)
    sig = torch.empty(B, device=device); rgb = torch.empty(B, 3, device=device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    out = {}

    def time_it(fn, iters=20):
        for _ in range(3):
            fn()
        evs = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b) for a, b in evs)
        return ts[len(ts) // 2] * 1e-3

    for name, xs, ds in (("random", x_rand, d), ("coherent", x_coh, d_coh)):
        t_f = time_it(lambda: field(xs, ds, out_sigmas=sig, out_rgbs=rgb))
        x01 = ((xs + 1) / 2).contiguous()
        feat = torch.empty(B, 32, dtype=torch.half, device=device)
        t_g = time_it(lambda: L.call("ntx_grid_encode_forward", L.ptr(x01), L.ptr(field.table), L.ptr(field.offsets), L.ptr(feat), B, 3, 2, 16, field.S,
                                     field.H, 0, None, 0, 1, L.F16, L.LAYOUT_BLC, L.stream()))
        out[name] = {"fused_field_msamples_per_s": B / t_f / 1e6, "fused_field_us": t_f * 1e6,
                     "fused_field_gbs": B * FIELD_BYTES_PER_SAMPLE / t_f / 1e9, "fused_field_frac_hbm": B * FIELD_BYTES_PER_SAMPLE / t_f / 1e9 / peaks["hbm_gbs"],
                     "fused_field_tflops": B * 36864 / t_f / 1e12,
                     "grid_encode_msamples_per_s": B / t_g / 1e6, "grid_encode_us": t_g * 1e6, "grid_encode_gbs": B * GRID_BYTES_PER_SAMPLE / t_g / 1e9,
                     "grid_encode_frac_hbm": B * GRID_BYTES_PER_SAMPLE / t_g / 1e9 / peaks["hbm_gbs"]}
    feat = torch.randn(B, 32, device=device).half()
    h = torch.empty(B, 16, dtype=torch.half, device=device)
    t_m = time_it(lambda: L.call("ntx_ffmlp_inference", L.ptr(feat), L.ptr(field.w_sigma), B, 32, 16, 64, 2, 0, 6, None, L.ptr(h), L.stream()))
    out["ffmlp_32_64_64_16"] = {"us": t_m * 1e6, "tflops": B * 14336 / t_m / 1e12, "frac_tensor_peak": B * 14336 / t_m / 1e12 / peaks["bf16_tflops"],
                                "io_gbs": B * 96 / t_m / 1e9, "io_frac_hbm": B * 96 / t_m / 1e9 / peaks["hbm_gbs"]}
    out["note"] = "2^20 samples, fp16 table 23.3 MiB (L2-resident), L2 flushed before every timed launch, median of 20"
    return out


if __name__ == "__main__":
    main()
