"""ctypes binding of the C-ABI library ``libnvsf_b200.so`` (include/nvsf_b200.h).

This is the whole "thin C-ABI torch-extension layer": tensors are passed as raw
device pointers plus the current CUDA stream handle; nothing torch-specific
crosses the boundary.  There is no fallback — if the library is missing or a
call fails the caller gets an exception.
"""
import ctypes
import contextlib
import functools
import threading
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# NVSF_B200_LIB: development override (A/B builds of the same sources); default = the in-tree library
LIB_PATH = os.environ.get("NVSF_B200_LIB") or os.path.join(_HERE, "libnvsf_b200.so")

_p = ctypes.c_void_p
_u32 = ctypes.c_uint32
_f32 = ctypes.c_float
_sz = ctypes.c_size_t
_int = ctypes.c_int

# name -> (restype, argtypes); mirrors include/nvsf_b200.h one to one.
PROTOTYPES = {
    "nvsf_abi_version": (_int, []),
    "nvsf_status_string": (ctypes.c_char_p, [_int]),
    "nvsf_near_far_from_aabb": (_int, [_p, _p, _p, _u32, _f32, _p, _p, _p]),
    "nvsf_sph_from_ray": (_int, [_p, _p, _f32, _u32, _p, _p]),
    "nvsf_morton3D": (_int, [_p, _u32, _p, _p]),
    "nvsf_morton3D_invert": (_int, [_p, _u32, _p, _p]),
    "nvsf_packbits": (_int, [_p, _u32, _f32, _p, _p]),
    "nvsf_march_rays_train_workspace_bytes": (_sz, [_u32]),
    "nvsf_march_rays_train": (
        _int,
        [_p, _p, _p, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _p, _p,
         _p, _sz, _p],
    ),
    "nvsf_march_rays_train_count": (
        _int,
        [_p, _p, _p, _f32, _f32, _u32, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _sz, _p],
    ),
    "nvsf_march_rays_train_write": (
        _int,
        [_p, _p, _p, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _p, _p,
         _u32, _p],
    ),
    "nvsf_march_rays_train_write_ws": (
        _int,
        [_p, _p, _p, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _p, _p,
         _u32, _p, _sz, _p],
    ),
    "nvsf_composite_rays_train_forward": (
        _int, [_p, _p, _p, _p, _u32, _u32, _f32, _p, _p, _p, _p]),
    "nvsf_composite_rays_train_backward": (
        _int, [_p, _p, _p, _p, _p, _p, _p, _p, _u32, _u32, _f32, _p, _p, _p]),
    "nvsf_march_rays": (
        _int,
        [_u32, _u32, _p, _p, _p, _p, _f32, _f32, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _p,
         _u32, _p],
    ),
    "nvsf_composite_rays": (_int, [_u32, _u32, _f32, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    # Part 2 (struct pointers are refined to typed pointers in field.py)
    "nvsf_field_workspace_bytes": (_sz, [_p]),
    "nvsf_field_pack_params": (_int, [_p, _p, _u32, _p, _sz, _p]),
    "nvsf_field_pack_time": (_int, [_p, _p, _p, _p, _sz, _p]),
    "nvsf_field_density_scratch_bytes": (_sz, [_u32]),
    "nvsf_field_density": (_int, [_p, _p, _p, _u32, _p, _p, _p, _p, _p, _sz, _p]),
    "nvsf_set_option": (_int, [ctypes.c_char_p, _int]),
    "nvsf_density_mode_get": (_int, []),
    "nvsf_get_option": (_int, [ctypes.c_char_p]),
    "nvsf_stage_timing_read": (_int, [_p, _p]),
    "nvsf_render_uniform_scratch_bytes": (_sz, [_u32, _u32]),
    "nvsf_render_uniform_density": (_int, [_p, _p, _p, _p, _p, _p, _p, _u32, _u32, _p, _sz, _p]),
    "nvsf_render_uniform_composite": (_int, [_p, _p, _u32, _p, _p, _p, _p, _u32, _u32, _f32, _p, _sz,
                                             _p, _p, _p, _p, _p, _p]),
    "nvsf_render_uniform": (_int, [_p, _p, _u32, _p, _p, _p, _p, _p, _u32, _u32, _f32, _p, _sz, _p,
                                   _p, _p, _p, _p, _p]),
    # Part 3 — training
    "nvsf_render_uniform_saved_bytes": (_sz, [_u32, _u32]),
    "nvsf_render_uniform_backward_scratch_bytes": (_sz, [_p, _u32, _u32]),
    "nvsf_render_uniform_debug_layout": (None, [_p, _u32, _u32, _p]),
    "nvsf_render_uniform_train_forward": (_int, [_p, _p, _u32, _p, _p, _p, _p, _p, _u32, _u32, _f32, _p,
                                                 _sz, _p, _p, _p, _p, _p, _p]),
    "nvsf_render_uniform_backward": (_int, [_p, _p, _p, _u32, _p, _p, _p, _p, _p, _u32, _u32, _f32, _p,
                                            _sz, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "nvsf_field_flow_scratch_bytes": (_sz, [_p, _u32]),
    "nvsf_field_flow_forward": (_int, [_p, _p, _p, _u32, _p, _p, _p, _sz, _p]),
    "nvsf_field_flow_backward": (_int, [_p, _p, _p, _p, _u32, _p, _p, _p, _p, _p, _sz, _p]),
    "nvsf_adam_step": (_int, [_p, _p, _p, _p, _sz, _f32, _f32, _f32, _f32, _u32, _f32, _p]),
    "nvsf_grad_found_inf": (_int, [_p, _sz, _p, _p]),
    "nvsf_adam_begin": (_int, [_p, _p, _f32, _f32, _p]),
    "nvsf_adam_step_guarded": (_int, [_p, _p, _p, _p, _sz, _f32, _f32, _f32, _f32, _p, _f32, _p]),
    "nvsf_ema_update": (_int, [_p, _p, _sz, _f32, _p]),
    "nvsf_field_color": (_int, [_p, _p, _u32, _p, _p, _u32, _u32, _p, _u32, _p, _u32, _p]),
    # Part 4 — ray generation, occupancy grid, alive-list compaction
    "nvsf_get_lidar_rays": (_int, [_p, _p, _u32, _u32, _u32, _f32, _f32, _f32, _p, _p, _p]),
    "nvsf_get_rays": (_int, [_p, _p, _u32, _u32, _u32, _f32, _f32, _f32, _f32, _p, _p, _p]),
    "nvsf_error_map_sample": (_int, [_p, _p, _p, _u32, _u32, _u32, _u32, _p, _p, _p]),
    "nvsf_error_map_update": (_int, [_p, _u32, _p, _u32, _p, _p]),
    "nvsf_grid_cell_points": (_int, [_u32, _u32, _f32, _p, _p, _p]),
    "nvsf_grid_cell_points_range": (_int, [_u32, _u32, _f32, _p, ctypes.c_uint64, ctypes.c_uint64, _p, _p]),
    "nvsf_grid_accumulate": (_int, [_p, _p, _u32, _f32, _u32, _p]),
    "nvsf_grid_update_workspace_bytes": (_sz, [_u32]),
    "nvsf_grid_update": (_int, [_p, _p, _u32, _f32, _f32, _p, _p, _p, _sz, _p]),
    "nvsf_compact_alive_workspace_bytes": (_sz, [_u32]),
    "nvsf_compact_alive": (_int, [_p, _u32, _p, _p, _p, _sz, _p]),
    # Part 5 — loss head
    "nvsf_loss_lidar": (_int, [_p, _p, _p, _u32, _p, _p, _p, _p, _p]),
    "nvsf_loss_elementwise": (_int, [_p, _p, _sz, _int, _f32, _f32, _p, _p, _p]),
    "nvsf_loss_los": (_int, [_p, _p, _p, _u32, _u32, _f32, _p, _p, _p, _sz, _p]),
    "nvsf_patch_grad_masks": (_int, [_p, _u32, _u32, _p, _u32, _u32, _u32, _f32, _f32, _p, _p, _p]),
    "nvsf_loss_patch": (_int, [_p, _p, _p, _p, _p, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _p]),
    "nvsf_chamfer_workspace_bytes": (_sz, [_u32, _u32, _u32]),
    "nvsf_chamfer_forward": (_int, [_p, _p, _u32, _u32, _u32, _p, _p, _p, _p, _p, _sz, _p]),
    "nvsf_chamfer_backward": (_int, [_p, _p, _u32, _u32, _u32, _p, _p, _p, _p, _p, _p, _p]),
    # Part 6 — evaluation
    "nvsf_chamfer_forward_counted": (_int, [_p, _p, _u32, _u32, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "nvsf_lidar_points_workspace_bytes": (_sz, [_u32, _u32]),
    "nvsf_lidar_points": (_int, [_p, _p, _f32, _p, _u32, _u32, _f32, _f32, _f32, _f32, _p, _p, _p, _sz, _p]),
    "nvsf_range_image_workspace_bytes": (_sz, [_u32, _u32, _u32]),
    "nvsf_range_image": (_int, [_p, _u32, _p, _u32, _u32, _p, _u32, _u32, _f32, _f32, _f32, _f32, _f32, _p, _p, _p,
                                _sz, _p]),
    "nvsf_eval_lidar_workspace_bytes": (_sz, [_u32, _u32]),
    "nvsf_eval_lidar": (_int, [_p, _p, _p, _u32, _u32, _f32, _f32, _f32, _f32, _f32, _f32, _p, _p, _sz, _p]),
    "nvsf_eval_camera_workspace_bytes": (_sz, [_u32, _u32]),
    "nvsf_eval_camera": (_int, [_p, _p, _u32, _u32, _p, _p, _sz, _p]),
    # Part 7 — mesh extraction
    "nvsf_marching_cubes_workspace_bytes": (_sz, [_u32, _u32, _u32]),
    "nvsf_marching_cubes_count": (_int, [_p, _u32, _u32, _u32, _f32, _p, _p, _sz, _p]),
    "nvsf_marching_cubes_write": (_int, [_p, _u32, _u32, _u32, _f32, _p, ctypes.c_uint64, _p, ctypes.c_uint64, _p,
                                         _sz, _p]),
}

_lib = None


class NvsfError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raise loudly if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA library has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`). "
            "nvsf_b200 has no CPU or PyTorch fallback."
        )
    handle = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(handle, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    got = handle.nvsf_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libnvsf_b200.so ABI {got} != python binding ABI {ABI_VERSION}; rebuild")
    _lib = handle
    return _lib


ABI_VERSION = 17


def check(status, what=""):
    if status != 0:
        msg = lib().nvsf_status_string(status).decode()
        raise NvsfError(f"{what}: {msg} (status {status})")


# ---- tuning options: process-wide in the C ABI, per model in this host mirror ----------------------------------
# nvsf_set_option writes process-wide switches that the launch code reads on the host at launch time.  The host
# mirror gives them per-model meaning and makes them safe with worker threads: every entry point of NeRFNetwork
# runs inside option_scope(model.options) — one re-entrant lock around "apply this model's overrides, enqueue the
# launches, restore" (the kernels themselves run asynchronously, outside the lock).
_OPTION_LOCK = threading.RLock()
_OPTION_LOCK_TIMEOUT_S = 120.0


def _acquire_option_lock():
    if not _OPTION_LOCK.acquire(timeout=_OPTION_LOCK_TIMEOUT_S):
        raise NvsfError(f"the option lock has been held by another thread for {_OPTION_LOCK_TIMEOUT_S:.0f} s "
                        "(is .backward() running inside a hand-opened option_scope? pass options=... to the model)")


@contextlib.contextmanager
def option_scope(overrides=None):
    """Hold the option lock; with `overrides` ({name: int}) set them for the duration and restore the previous
    values afterwards.  Unknown names / rejected values raise NvsfError before anything is launched."""
    # (a bounded wait: a thread that opens a scope by hand and calls loss.backward() inside it would otherwise wait
    #  forever for the autograd thread, which needs the same lock — give the MODEL its options instead)
    _acquire_option_lock()
    try:
        if not overrides:
            yield
            return
        L = lib()
        saved = []
        try:
            for name, value in overrides.items():
                key = name.encode()
                old = L.nvsf_get_option(key)
                check(L.nvsf_set_option(key, int(value)), f"set_option({name}={value})")
                saved.append((key, old))
            yield
        finally:
            for key, old in reversed(saved):
                L.nvsf_set_option(key, old)
    finally:
        _OPTION_LOCK.release()


def with_options(fn):
    """Method decorator: run under option_scope(self.options) (see above)."""

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with option_scope(getattr(self, "options", None)):
            return fn(self, *args, **kwargs)

    return wrapper


def ptr(t):
    """Raw device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr() or None


def stream_ptr():
    import torch

    return torch.cuda.current_stream().cuda_stream or None


def device_guard(fn):
    """Run `fn` with the CUDA device of its first CUDA tensor (or of the first nn.Module with CUDA
    parameters) current, as torch's own extensions do through their device guard: the kernels behind
    the C ABI launch on the current device and on its current stream (`stream_ptr`)."""
    import torch

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        for a in args:
            if isinstance(a, torch.Tensor):
                if a.is_cuda:
                    dev = a.device
                    break
            elif isinstance(a, torch.nn.Module):
                p = next(a.parameters(), None)
                if p is not None and p.is_cuda:
                    dev = p.device
                    break
        # the option lock: a launch never observes another thread's model-scoped overrides half applied
        _acquire_option_lock()
        try:
            if dev is None or dev.index == torch.cuda.current_device():
                return fn(*args, **kwargs)
            with torch.cuda.device(dev):
                return fn(*args, **kwargs)
        finally:
            _OPTION_LOCK.release()

    return wrapper
