"""ctypes binding of libntx.so (the C ABI declared in include/ntx.h).

There is deliberately no CPU fallback: if the library is missing or a call fails, a RuntimeError is raised —
the same exception type the reference's TORCH_CHECK / std::runtime_error surface as in Python.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NTX_LIB_PATH") or os.path.join(_HERE, "lib", "libntx.so")   # NTX_LIB_PATH: development (tools/tune.py variants)
_lib = None

F32, F16, F64 = 0, 1, 2
LAYOUT_LBC, LAYOUT_BLC = 0, 1
_DTYPE_ID = {torch.float32: F32, torch.float16: F16, torch.float64: F64}

_u32, _f32, _int, _vp, _sz = C.c_uint32, C.c_float, C.c_int, C.c_void_p, C.c_size_t
_SIGS = {
    "ntx_grid_encode_forward": [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _f32, _u32, _int, _vp, _u32, _int, _int, _int, _vp],
    "ntx_grid_encode_backward": [_vp, _vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _f32, _u32, _int, _vp, _vp, _u32, _int, _int, _int, _vp],
    "ntx_grid_level_scales": [_f32, _u32, _u32, _vp, _vp],
    "ntx_grid_debug_indices": [_vp, _vp, _u32, _u32, _u32, _f32, _u32, _u32, _int, _vp, _vp],
    "ntx_ffmlp_forward": [_vp, _vp, _u32, _u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp],
    "ntx_ffmlp_inference": [_vp, _vp, _u32, _u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp],
    "ntx_ffmlp_backward": [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _u32, _u32, _u32, _int, _vp, _vp, _vp, _vp, _vp],
    "ntx_allocate_splitk": [_sz],
    "ntx_free_splitk": [],
    "ntx_sh_encode_forward": [_vp, _vp, _u32, _u32, _u32, _int, _vp, _vp],
    "ntx_sh_encode_backward": [_vp, _vp, _u32, _u32, _u32, _vp, _vp, _vp],
    "ntx_near_far_from_aabb": [_vp, _vp, _vp, _u32, _f32, _vp, _vp, _vp],
    "ntx_polar_from_ray": [_vp, _vp, _f32, _u32, _vp, _vp],
    "ntx_morton3D": [_vp, _u32, _vp, _vp],
    "ntx_morton3D_invert": [_vp, _u32, _vp, _vp],
    "ntx_packbits": [_vp, _u32, _f32, _vp, _vp],
    "ntx_march_rays_train": [_vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _vp, _vp],
    "ntx_composite_rays_train_forward": [_vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp],
    "ntx_composite_rays_train_backward": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp],
    "ntx_march_rays": [_u32, _u32, _vp, _vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _int, _u32, _vp, _vp],
    "ntx_build_occupancy_mip": [_vp, _u32, _u32, _vp, _vp],
    "ntx_composite_rays": [_u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "ntx_compact_rays": [_u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "ntx_ngp_field_forward": [_vp, _vp, _vp, _u32, _f32, _vp, _vp, _u32, _f32, _u32, _int, _vp, _vp, _f32, _vp, _vp, _vp],
    "ntx_render_rays": [_vp, _vp, _u32, _vp, _f32, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _u32, _f32, _u32, _int, _vp, _vp, _f32,
                        _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "ntx_unshard_frame": [_vp, _u32, _u32, _u32, _u32, _f32, _vp, _vp, _vp, _vp],
    "ntx_unshard_frame_peers": [_vp, _sz, _u32, _u32, _u32, _u32, _f32, _vp, _vp, _vp, _vp],
    "ntx_mesh_create": [_vp, _u32, _vp, _u32, _vp],
    "ntx_mesh_destroy": [_vp],
    "ntx_mesh_info": [_vp, _vp],
    "ntx_mesh_trace": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _vp],
    "ntx_mesh_knn": [_vp, _vp, _u32, _u32, _f32, _vp, _vp, _vp],
    "ntx_mesh_project": [_vp, _vp, _vp, _u32, _u32, _f32, _f32, _vp, _vp, _vp, _vp, _vp],
    "ntx_texture_field_density": [_vp, _vp, _vp, _u32, _u32, _f32, _f32, _f32, _f32, _vp, _vp, _u32, _f32, _u32, _int, _vp, _vp, _vp, _vp],
    "ntx_update_density_grid": [_vp, _vp, _u32, _u32, _f32, _f32, _f32, _f32, _vp, _vp, _u32, _f32, _u32, _int, _vp, _vp, _u32, _vp, _int, _vp, _vp, _vp],
}
_SIZE_FNS = {
    "ntx_update_density_grid_workspace_bytes": [_u32, _u32],
    "ntx_march_rays_train_workspace_bytes": [_u32],
    "ntx_compact_rays_workspace_bytes": [_u32],
    "ntx_occupancy_mip_bytes": [_u32, _u32],
    "ntx_render_rays_workspace_bytes": [_u32, _u32],
    "ntx_ffmlp_backward_workspace_bytes": [_u32, _u32, _u32, _u32],
}


def lib():
    """Load libntx.so (building is the job of __graft_entry__.build() / `python -m nerf_texture_b200.build`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libntx.so not found at %s — build it with `python -m nerf_texture_b200.build` (there is no CPU fallback)" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        l.ntx_last_error.restype = C.c_char_p
        for name, sig in _SIGS.items():
            if hasattr(l, name):
                fn = getattr(l, name)
                fn.argtypes = sig
                fn.restype = C.c_int
        for name, sig in _SIZE_FNS.items():
            if hasattr(l, name):
                fn = getattr(l, name)
                fn.argtypes = sig
                fn.restype = C.c_size_t
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError(lib().ntx_last_error().decode() or "libntx error %d" % rc)


launches = 0  # number of libntx kernel-launching calls made by this process (bench.py reports the delta as gpu_launches)
_NO_LAUNCH = {"ntx_allocate_splitk", "ntx_free_splitk", "ntx_mesh_create", "ntx_mesh_destroy", "ntx_mesh_info"}


def call(name, *args):
    global launches
    check(getattr(lib(), name)(*args))
    if name not in _NO_LAUNCH:
        launches += 1


def ptr(t, dtype=None):
    """device pointer of a CUDA tensor (None -> NULL); the reference's CHECK_CUDA / CHECK_CONTIGUOUS / CHECK_IS_INT /
    CHECK_IS_FLOATING live here: a wrong dtype or a tensor on another GPU raises instead of being reinterpreted
    (the reference raises through data_ptr<T>() in that case)"""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("tensor must be a CUDA tensor")
    if not t.is_contiguous():
        raise RuntimeError("tensor must be a contiguous tensor")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("tensor must be a %s tensor (got %s)" % (str(dtype).replace("torch.", ""), str(t.dtype).replace("torch.", "")))
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError("tensor is on cuda:%d but the current device is cuda:%d" % (t.device.index, torch.cuda.current_device()))
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def dtype_id(dt):
    if dt not in _DTYPE_ID:
        raise RuntimeError("tensor must be a floating tensor")
    return _DTYPE_ID[dt]


_workspaces = {}


def workspace(kind, nbytes, device):
    """Zero-initialised, self-cleaning scan workspace, one per (kind, device, stream) and grown on demand."""
    key = (kind, device.index, stream())
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(int(nbytes), 4096), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def bind_host_thread_to_gpu(device_index):
    """Pin the calling thread (and what it allocates next: pinned staging buffers, the frame mailbox) to the CPUs of the NUMA node the
    GPU hangs off (NVML's ideal CPU affinity).  On a two-socket B200 box a rank whose pinned buffers live on the far socket pays for it
    in every host<->device copy and every mailbox read; returns the previous affinity (for os.sched_setaffinity) or None if NVML is
    not available.  Best effort: never raises."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        prev = os.sched_getaffinity(0)
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(int(device_index)))
        return prev
    except Exception:
        return None
