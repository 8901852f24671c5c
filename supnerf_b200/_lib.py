"""ctypes binding of libsupnerf_b200.so (the C ABI declared in include/supnerf_b200.h).

There is no fallback: if the library is missing, or a call fails, this raises."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsupnerf_b200.so")

c_f = ctypes.c_void_p  # device float*
c_i64, c_i32, c_flt, c_sz = ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_size_t


class SnbArch(ctypes.Structure):
    _fields_ = [("arch", c_i32), ("shape_blocks", c_i32), ("texture_blocks", c_i32), ("W", c_i32),
                ("latent_dim", c_i32), ("num_xyz_freq", c_i32), ("num_dir_freq", c_i32)]


class SnbRenderDesc(ctypes.Structure):
    _fields_ = [("n_rays", c_i64), ("n_samples", c_i32), ("precision", c_i32), ("flags", c_i32), ("half_diag", c_flt),
                ("aabb_half", c_flt * 3), ("mode", c_i32), ("obj_diag", c_flt), ("shapenet_swap", c_i32)]


class SnbBatchDesc(ctypes.Structure):
    _fields_ = [("n_objs", c_i32), ("n_samples", c_i32), ("rays_per_obj", c_i64), ("flags", c_i32), ("reserved", c_i32)]


class SnbShellBatchDesc(ctypes.Structure):
    _fields_ = [("n_objs", c_i32), ("n_samples", c_i32), ("rays_per_obj", c_i64), ("precision", c_i32), ("flags", c_i32),
                ("shapenet_swap", c_i32), ("reserved", c_i32)]


# name -> (restype, argtypes); mirrors include/supnerf_b200.h one to one
SIGNATURES = {
    "snb_abi_version": (c_i32, []),
    "snb_last_error": (ctypes.c_char_p, []),
    "snb_launch_count": (ctypes.c_uint64, []),
    "snb_device_info": (c_i32, [ctypes.POINTER(c_i32)] * 3),
    "snb_composite_fwd": (c_i32, [c_f, c_f, c_f, c_i64, c_i64, c_i32, c_i32, c_f, c_f, c_f, c_f]),
    "snb_composite_bwd": (c_i32, [c_f, c_f, c_f, c_i64, c_i64, c_i32, c_i32, c_f, c_f, c_f, c_f, c_f, c_f, c_f]),
    "snb_get_rays_fwd": (c_i32, [c_f, c_f, c_i64, c_f, c_f, c_f, c_f, c_f]),
    "snb_get_rays_bwd": (c_i32, [c_f, c_f, c_i64, c_f, c_f, c_f, c_f, c_f, c_f]),
    "snb_ray_box_fwd": (c_i32, [c_f, c_f, c_f, c_f, c_i64, c_f, c_f, c_f, c_f]),
    "snb_ray_box_bwd": (c_i32, [c_f, c_f, c_f, c_f, c_i64, c_f, c_f, c_f, c_f, c_f, c_f, c_f]),
    "snb_sample_box_fwd": (c_i32, [c_f, c_f, c_f, c_f, c_i64, c_i32, c_flt, ctypes.POINTER(c_flt), c_f, c_f, c_f, c_f, c_f]),
    "snb_sample_box_bwd": (c_i32, [c_f, c_f, c_f, c_f, c_i64, c_i32, c_flt, ctypes.POINTER(c_flt), c_f, c_f, c_f, c_f, c_f, c_i32, c_f]),
    "snb_stratified_z_fwd": (c_i32, [c_f, c_i32, c_f, c_f, c_i64, c_i32, c_f, c_f]),
    "snb_stratified_z_bwd": (c_i32, [c_f, c_f, c_i64, c_i32, c_f, c_f, c_f, c_f]),
    "snb_sample_shell_fwd": (c_i32, [c_f, c_f, c_f, c_i64, c_i32, c_flt, c_i32, c_f, c_f, c_f]),
    "snb_sample_shell_bwd": (c_i32, [c_f, c_i64, c_i32, c_flt, c_i32, c_f, c_f, c_f, c_f, c_f]),
    "snb_jitter_fill": (c_i32, [ctypes.c_uint64, c_f, c_i64, c_i32, c_f, c_f]),
    "snb_create": (c_i32, [ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(SnbArch)]),
    "snb_destroy": (c_i32, [ctypes.c_void_p]),
    "snb_num_weight_tensors": (c_i32, [ctypes.c_void_p]),
    "snb_layer_shape": (c_i32, [ctypes.c_void_p, c_i32, ctypes.POINTER(c_i32), ctypes.POINTER(c_i32)]),
    "snb_set_weights": (c_i32, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), c_i32]),
    "snb_packed_bytes": (c_sz, [ctypes.c_void_p]),
    "snb_tc_set_debug": (c_i32, [ctypes.c_void_p, c_f]),
    "snb_tc_set_trace": (c_i32, [ctypes.c_void_p, c_f]),
    "snb_tc_set_cg2": (c_i32, [ctypes.c_void_p, c_i32]),
    "snb_kernel_timing_enable": (c_i32, [ctypes.c_void_p, c_i32]),
    "snb_kernel_timing_read": (c_i32, [ctypes.c_void_p, c_i32, ctypes.POINTER(c_flt), c_i32]),
    "snb_pack_weights": (c_i32, [ctypes.c_void_p, c_f, c_f]),
    "snb_mlp_workspace_bytes": (c_sz, [ctypes.c_void_p, c_i64, c_i64, c_i32]),
    "snb_mlp_bwd_scratch_bytes": (c_sz, [ctypes.c_void_p, c_i64, c_i64, c_i32]),
    "snb_mlp_fwd": (c_i32, [ctypes.c_void_p, c_i32, c_f, c_f, c_i64, c_i64, c_f, c_f, c_f, c_f, c_f, c_f]),
    "snb_mlp_bwd": (c_i32, [ctypes.c_void_p, c_i32, c_f, c_f, c_i64, c_i64, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_f,
                            c_f, c_f, ctypes.POINTER(ctypes.c_void_p), c_f]),
    "snb_refine_loss_scratch_bytes": (c_sz, []),
    "snb_refine_loss_fwd": (c_i32, [c_f, c_f, c_f, c_f, c_i64, c_flt, c_f, c_f, c_f, c_f]),
    "snb_refine_loss_bwd": (c_i32, [c_f, c_f, c_f, c_f, c_i64, c_flt, c_f, c_f, c_f, c_f, c_f]),
    "snb_merge_sort_samples": (c_i32, [c_f, c_f, c_f, c_i64, c_i32, c_f, c_f, c_f, c_f, c_f]),
    "snb_render_workspace_bytes": (c_sz, [ctypes.c_void_p, ctypes.POINTER(SnbRenderDesc)]),
    "snb_render_bwd_scratch_bytes": (c_sz, [ctypes.c_void_p, ctypes.POINTER(SnbRenderDesc)]),
    "snb_render_fwd": (c_i32, [ctypes.c_void_p, ctypes.POINTER(SnbRenderDesc)] + [c_f] * 14),
    "snb_render_bwd": (c_i32, [ctypes.c_void_p, ctypes.POINTER(SnbRenderDesc)] + [c_f] * 16 + [ctypes.POINTER(ctypes.c_void_p), c_f]),
    "snb_allreduce_grads": (c_i32, [ctypes.c_void_p, ctypes.c_void_p, c_f, c_sz, c_f]),
    "snb_render_batch_workspace_bytes": (c_sz, [ctypes.c_void_p, ctypes.POINTER(SnbBatchDesc)]),
    "snb_render_batch_scratch_bytes": (c_sz, [ctypes.c_void_p, ctypes.POINTER(SnbBatchDesc)]),
    "snb_render_batch_fwd": (c_i32, [ctypes.c_void_p, ctypes.POINTER(SnbBatchDesc)] + [c_f] * 15),
    "snb_render_batch_bwd": (c_i32, [ctypes.c_void_p, ctypes.POINTER(SnbBatchDesc)] + [c_f] * 18),
    "snb_prepare_samples_batch": (c_i32, [c_f, c_f, c_f, c_f, c_f, c_f, c_f, c_i32, c_i64, c_i32, c_i32, c_f, c_f, c_f]),
    "snb_refine_loss_batch_scratch_bytes": (c_sz, [c_i32]),
    "snb_refine_loss_batch_fwd": (c_i32, [c_f, c_f, c_f, c_f, c_i32, c_i64, c_flt, c_f, c_f, c_f]),
    "snb_refine_loss_batch_bwd": (c_i32, [c_f, c_f, c_f, c_f, c_i32, c_i64, c_flt, c_f, c_f, c_f, c_f, c_f]),
    "snb_refine_pose_batch_bwd": (c_i32, [c_f, c_f, c_i32, c_i32, c_f, c_f, c_f, c_f]),
    "snb_refine_pose_slots_fwd": (c_i32, [c_f, c_f, c_i32, c_i32, c_f, c_i32, c_f, c_f, c_f, c_i32, c_f, c_f, c_f, c_f, c_f, c_f]),
    "snb_adamw_step_rows": (c_i32, [c_i32, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                    ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(c_i32), ctypes.POINTER(c_flt), c_flt, c_flt, c_flt, c_flt,
                                    c_i32, c_f, c_f, c_f, c_f, c_i32, c_f, c_i32, c_f]),
    "snb_render_shell_batch_workspace_bytes": (c_sz, [ctypes.c_void_p, ctypes.POINTER(SnbShellBatchDesc)]),
    "snb_render_shell_batch_scratch_bytes": (c_sz, [ctypes.c_void_p, ctypes.POINTER(SnbShellBatchDesc)]),
    "snb_render_shell_batch_fwd": (c_i32, [ctypes.c_void_p, ctypes.POINTER(SnbShellBatchDesc)] + [c_f] * 13),
    "snb_render_shell_batch_bwd": (c_i32, [ctypes.c_void_p, ctypes.POINTER(SnbShellBatchDesc)] + [c_f] * 17),
}

_lib = None


def load():
    """Load the shared library (once).  Raises if it has not been built — there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m supnerf_b200.build` (or __graft_entry__.build()). "
            "supnerf_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.snb_abi_version() != 2:
        raise ImportError("libsupnerf_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


class SnbError(RuntimeError):
    pass


def check(rc, what):
    if rc != 0:
        raise SnbError(f"{what} failed (rc={rc}): {load().snb_last_error().decode(errors='replace')}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  Tensors must be CUDA, fp32/uint8, contiguous."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    """cudaStream_t of torch's current stream on the current device (the raw accessor: torch.cuda.current_stream() builds a
    Stream object per call, ~10x the cost, and every C-ABI call needs this)."""
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NO_GUARD = _NoGuard()


def on_device(dev):
    """`with on_device(t.device):` == `with torch.cuda.device(t.device):`, but free when that device is already current."""
    if dev.index is None or torch._C._cuda_getDevice() == dev.index:
        return _NO_GUARD
    return torch.cuda.device(dev)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise SnbError("supnerf_b200 kernels need CUDA tensors; there is no CPU fallback")


def f32c(t):
    """contiguous fp32 view/copy on the same device"""
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()
