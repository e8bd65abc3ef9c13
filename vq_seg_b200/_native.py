"""ctypes binding of libvqseg.so (C ABI declared in include/vqseg.h).

There is NO CPU fallback: if the shared library is missing or the device is not a B200 the
calls raise.  Build with `python -m vq_seg_b200.build` (or `__graft_entry__.build()`).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvqseg.so")
DEV_LIB_PATH = os.path.join(_HERE, "libvqseg_dev.so")      # developer build (-DVQSEG_DEV): pipeline trace hooks, never shipped
_lib = None

i64, f32, vp, sz, ci = ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int

# name -> (restype, argtypes); mirrors include/vqseg.h one to one
SIGNATURES = {
    "vqseg_version": (ci, []),
    "vqseg_error_string": (ctypes.c_char_p, [ci]),
    "vqseg_codebook_blob_bytes": (sz, [i64, i64]),
    "vqseg_codebook_prepare_f32": (ci, [vp, i64, i64, vp, sz, vp]),
    "vqseg_codebook_prepare_ip_f32": (ci, [vp, i64, i64, vp, sz, vp]),
    "vqseg_samples_blob_bytes": (sz, [i64, i64]),
    "vqseg_samples_prepare_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, sz, vp]),
    "vqseg_assign_prepared_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, vp, i64, vp, vp, vp, ci, vp, sz, vp, vp]),
    "vqseg_assign_workspace_bytes": (sz, [i64, i64, i64, ci]),
    "vqseg_assign_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, vp, vp, vp, vp, i64, ci, ci, vp, sz, vp, vp]),
    "vqseg_unpack_keys": (ci, [vp, i64, vp, vp, vp, i64, vp]),
    "vqseg_gather_workspace_bytes": (sz, [i64, i64]),
    "vqseg_gather_ste_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, vp, vp, i64, i64, i64, vp, ci, vp, sz, vp]),
    "vqseg_forward_workspace_bytes": (sz, [i64, i64, i64]),
    "vqseg_vq_forward_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, vp, vp, vp, vp, vp, i64, i64, i64, vp,
                                  ci, ci, ci, vp, sz, vp, vp]),
    "vqseg_ste_bwd_f32": (ci, [vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64, vp, f32,
                               vp, i64, i64, i64, i64, i64, i64, vp]),
    "vqseg_rotate_bwd_f32": (ci, [vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64, vp, f32,
                                  vp, i64, i64, i64, i64, i64, i64, vp]),
    "vqseg_gather_bwd_codebook_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, vp, i64, vp]),
    "vqseg_code_stats_workspace_bytes": (sz, [i64, i64, i64, ci]),
    "vqseg_code_stats_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, vp, vp, ci, vp, sz, vp]),
    "vqseg_kmeans_finalize_f32": (ci, [vp, vp, vp, i64, i64, ci, vp]),
    "vqseg_code_usage": (ci, [vp, i64, vp, vp]),
    "vqseg_gather_rows_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, vp, vp]),
    "vqseg_l2norm_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, i64, i64, vp]),
    "vqseg_ema_update_f32": (ci, [vp, vp, vp, vp, vp, i64, i64, f32, f32, vp, vp]),
    "vqseg_ema_expire_workspace_bytes": (sz, [i64]),
    "vqseg_ema_update_expire_f32": (ci, [vp, vp, vp, vp, vp, i64, i64, f32, f32, f32, f32, vp, vp, vp, sz, vp]),
    "vqseg_dist_map_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, ci, vp, i64, i64, i64, vp, vp, vp, vp]),
    "vqseg_dist_map_bwd_f32": (ci, [vp, vp, i64, i64, i64, vp, i64, i64, i64, i64, i64, i64, vp, i64,
                                    vp, i64, i64, i64, vp, vp, vp]),
    "vqseg_sim_map_bwd_f32": (ci, [vp, i64, i64, i64, vp, i64, i64, i64, i64, i64, i64, vp, i64, vp, i64, i64, i64, vp, vp]),
    "vqseg_seghead_map_f32": (ci, [vp, i64, i64, i64, i64, i64, i64, vp, i64, ci, vp, i64, i64, i64, vp, vp, vp, ci, vp]),
    "vqseg_seghead_map_bwd_workspace_bytes": (sz, [i64, i64, i64, ci]),
    "vqseg_seghead_map_bwd_f32": (ci, [vp, vp, i64, i64, i64, vp, i64, i64, i64, i64, i64, i64, vp, i64, ci, vp,
                                       vp, i64, i64, i64, vp, ci, vp, sz, vp]),
}


class NativeLibraryError(RuntimeError):
    pass


def lib():
    """Loads libvqseg.so once; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                f"{LIB_PATH} not found: build it with `python -m vq_seg_b200.build`. "
                "vq_seg_b200 has no CPU / PyTorch fallback for its kernels.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError if the .so does not export it
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def use_dev_library():
    """scripts/gpu_dev.py only: bind the developer build (same ABI + vqseg_debug_set_trace) instead of the product .so."""
    global _lib
    handle = ctypes.CDLL(DEV_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)
        fn.restype, fn.argtypes = res, args
    handle.vqseg_debug_set_trace.restype, handle.vqseg_debug_set_trace.argtypes = None, [vp]
    _lib = handle
    return handle


class ProfileEvents:
    """Four caller-owned CUDA events handed to vqseg_assign_f32 / vqseg_vq_forward_f32 (`prof_events`): the call
    records [0],[1] around the tensor-core filter kernel and [2],[3] around the rescoring kernel."""

    def __init__(self):
        import torch
        self.events = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        for e in self.events:
            e.record()                      # torch creates the cudaEvent_t lazily, on the first record
        torch.cuda.synchronize()
        self.array = (vp * 4)(*[e.cuda_event for e in self.events])

    def _ms(self, a, b):
        try:                                # the caller has synchronised the stream / device
            return self.events[a].elapsed_time(self.events[b])
        except RuntimeError:
            return -1.0

    def filter_ms(self):
        return self._ms(0, 1)

    def rescore_ms(self):
        return self._ms(2, 3)


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().vqseg_error_string(rc).decode()
        raise RuntimeError(f"libvqseg {what} failed ({rc}): {msg}")
