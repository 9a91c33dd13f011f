"""Builds nerf_texture_b200/lib/libntx.so — the C-ABI CUDA library — with nvcc for sm_100a, in-tree.

    python -m nerf_texture_b200.build [--force] [--verbose]

Each .cu is compiled to an object (in parallel) and linked into one shared library with a static cudart, so the
.so only needs the CUDA driver on the GPU box.  No torch headers are involved: the kernels take raw pointers.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
# development variants: NTX_BUILD_TAG=probe NTX_NVCC_EXTRA=-DNTX_DEV_PROBES builds lib/libntx_probe.so next to the product library
# (select it at run time with NTX_LIB_PATH); the product build has no tag
_TAG = os.environ.get("NTX_BUILD_TAG", "")
OBJDIR = os.path.join(LIBDIR, "obj" + ("_" + _TAG if _TAG else ""))
LIB = os.path.join(LIBDIR, "libntx" + ("_" + _TAG if _TAG else "") + ".so")
# longest compile first (mlp.cu: ~55 s of ~100 s in all), so that a build with fewer jobs than sources is not left waiting on it at the end
SOURCES = ["mlp.cu", "grid.cu", "mlp_bwd.cu", "mesh.cu", "texture_field.cu", "raymarch.cu", "field.cu", "sh.cu", "api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr", "-Xptxas", "-v",
] + os.environ.get("NTX_NVCC_EXTRA", "").split()   # development only, e.g. -DNTX_DEV_PROBES (tools/field_probe.py)


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _deps(src):
    deps = [os.path.join(CSRC, src), os.path.join(HERE, "..", "include", "ntx.h")]
    deps += [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))]
    return deps


def _stamp(src):
    h = hashlib.sha1(" ".join(NVCC_FLAGS).encode())
    for d in sorted(_deps(src)):
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _compile(src, force, verbose):
    obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
    stamp_file = obj + ".stamp"
    stamp = _stamp(src)
    if not force and os.path.exists(obj) and os.path.exists(stamp_file) and open(stamp_file).read() == stamp:
        return obj, False, ""
    cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout[-6000:], r.stderr[-12000:]))
    with open(stamp_file, "w") as f:
        f.write(stamp)
    with open(obj + ".ptxas.log", "w") as f:
        f.write(r.stderr)
    return obj, True, r.stderr


def _mem_available_bytes():
    """memory this process can still use: MemAvailable, or less under a cgroup (v2) memory limit; None if unknown"""
    avail = None
    try:
        with open("/proc/meminfo") as f:
            avail = next(int(l.split()[1]) * 1024 for l in f if l.startswith("MemAvailable:"))
    except (OSError, StopIteration, ValueError):
        pass
    try:
        with open("/sys/fs/cgroup/memory.max") as f:
            limit = f.read().strip()
        if limit != "max":
            with open("/sys/fs/cgroup/memory.current") as f:
                free = int(limit) - int(f.read().strip())
            avail = free if avail is None else min(avail, free)
    except (OSError, ValueError):
        pass
    return avail


def _jobs(n):
    """parallel nvcc jobs: no more than the CPUs this process may run on (os.cpu_count() counts the host's in a container) and one per
    GB of available memory (cicc + ptxas of mlp.cu peak at ~0.6 GB, the other sources at ~0.25 GB)"""
    try:
        cpus = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        cpus = os.cpu_count() or 4
    mem = _mem_available_bytes()
    by_mem = max(1, mem // (1 << 30)) if mem is not None else cpus
    return max(1, min(n, cpus, by_mem))


def build(force=False, verbose=False):
    os.makedirs(OBJDIR, exist_ok=True)
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    with ThreadPoolExecutor(max_workers=_jobs(len(srcs))) as ex:
        results = list(ex.map(lambda s: _compile(s, force, verbose), srcs))
    objs = [r[0] for r in results]
    rebuilt = any(r[1] for r in results)
    if verbose:
        for s, r in zip(srcs, results):
            if r[1]:
                print("== %s ==\n%s" % (s, r[2]))
    if rebuilt or not os.path.exists(LIB):
        cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-cudart", "static", "-Xcompiler", "-fPIC"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv or "-v" in sys.argv))
